"""Read sets planned against the slot index's own geometry, so that its probe walks reach their edges on purpose.

TEST INFRASTRUCTURE.  Every stage reaches the prefix/suffix table through an open-addressing walk over 4-slot sectors that
starts in the key's home sector, moves on while a sector is full and wraps from the last sector of the index (or of the
key's shard) to its first.  A random key homes in the last sector with probability 1 / nsec, so the ordinary data sets wrap
and build long chains only by chance.  The sets here fix the number of unique reads U first, which fixes the index size
(table_shard_slots in csrc/table.cu, restated below), and then choose keys by rejection sampling so that they home where a
chain has to form:

  wrap_end      the last 8 sectors of the single table overfilled: the chain runs past nsec - 1 and on from sector 0
  long_run      16 or more consecutive full sectors in the middle of the index: one read probes a long walk and short ones
  bucket_seam   a chain across the boundary between two slot ranges of the bucketed build (a bucket = top 8 hash bits)
  shard_ends2/3 chains that wrap at the end of shard 0 and of shard 1 of a 2- / 3-shard table

Hashes, home sectors, owners and tags come from tests/table_ref.py, which restates core.cuh.

The crafted keys sit in a genome: block j of D bases is the crafted h-mer (or its reverse complement) and a random spacer.
The read of block j starts at the block (forward) or ends at its h-mer (a reverse-strand read, given reverse complemented),
and two spacer bases are fixed to A so that every crafted read is stored in the orientation planned: its first h bases are
then the key of the type planned (0 / 2 as given, 1 / 3 through their reverse complement).  A read spans the next block's
h-mer too, and a second read starts 7 bases into every block, so the crafted keys are also interior windows of the search.
A masked key (110 reads) and a run key (40 reads) share their first h bases with distinct remainders and home at the end of
the crowded chain with the largest hashes of their sector, so that the reference build (keys in hash order) puts them in
the part of the chain that was pushed furthest (past the wrap where there is one).  Random reads fill the set up to U.
"""
from __future__ import annotations

import functools

import numpy as np

import table_ref

SETS = ["wrap_end", "long_run", "bucket_seam", "shard_ends2", "shard_ends3"]
KS = [32, 45, 70]
U_PLAN = 3000
MASKED_READS, RUN_READS = 110, 40
BUCKET = 128                         # bucket_seam: the chain crosses from bucket 127 into bucket 128
LONG_RUN_SECTORS, LONG_WALK = 16, 10
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_u = np.uint64

# (block length D, read length L) per h: the last base of a forward read and the first base of a reverse-strand read fall in
# the spacer of a block ((L - 1) % D and (h - L) % D are both >= h), and a read spans the next block's h-mer (D + h <= L)
GEOMETRY = {32: (50, 100), 45: (60, 120), 64: (80, 150)}


def table_sectors(U: int, world: int = 1) -> int:
    """sectors of one shard of the slot index (csrc/table.cu table_shard_slots)"""
    n = 4 * U
    nsec = (n + n // 2 + 3) // 4
    if world > 1:
        nsec = nsec // world + nsec // (10 * world) + 1
    return max(nsec, 256)


def world_of(name: str) -> int:
    return int(name[-1]) if name.startswith("shard_ends") else 1


def _key_words(codes: np.ndarray, h: int):
    """(v0, v1) of h-mers given as rows of 2-bit codes (table_ref.Keys' fold)"""
    w = codes.astype(np.uint64)
    v0 = np.zeros(len(codes), np.uint64)
    v1 = np.zeros(len(codes), np.uint64)
    split = max(h - 32, 0)
    for t in range(split):
        v0 = (v0 << _u(2)) | w[:, t]
    for t in range(split, h):
        v1 = (v1 << _u(2)) | w[:, t]
    return v0, v1


def _hash(codes: np.ndarray, h: int) -> np.ndarray:
    return table_ref.hash_key(*_key_words(codes, h))


def _rc(codes: np.ndarray) -> np.ndarray:
    return (3 - codes)[..., ::-1]


class _Sampler:
    """h-mers drawn in batches of random candidates; a draw takes the first unused candidate that meets its target"""

    def __init__(self, rng, h, nsec, world):
        self.rng, self.h, self.nsec, self.world = rng, h, nsec, world
        self.pools = {}

    def _pool(self, first, target_rc):
        if (first, target_rc) not in self.pools:
            c = self.rng.integers(0, 4, size=(400_000, self.h), dtype=np.uint8)
            c[:, 0] = first
            hsh = _hash(_rc(c) if target_rc else c, self.h)
            with np.errstate(over="ignore"):      # an eighth of a sector further is the next sector (or past 2^64)
                up = hsh + _u(1 << 61) // _u(self.nsec)
            sec = table_ref.home_sector(hsh, self.nsec).astype(np.int64)
            top = (up < hsh) | (table_ref.home_sector(up, self.nsec).astype(np.int64) > sec)
            self.pools[first, target_rc] = [c, hsh, sec, top, table_ref.key_owner(hsh, self.world), np.zeros(len(c), bool)]
        return self.pools[first, target_rc]

    def draw(self, first: int, target_rc: bool, lo: int, hi: int, owner: int = 0, top: bool = False):
        """an h-mer starting with base `first` whose key (its reverse complement when target_rc) homes in [lo, hi) of the
        shard `owner`; top: in the top eighth of its home sector's hash range"""
        c, hsh, sec, is_top, own, used = self._pool(first, target_rc)
        ok = (sec >= lo) & (sec < hi) & (own == owner) & ~used
        if top:
            ok &= is_top
        at = np.flatnonzero(ok)
        assert len(at), "no h-mer found for the target"
        used[at[0]] = True
        return c[at[0]]


class Plan:
    """A planned set: reads (bytes, as given to the pipeline), k, h, U, world, nsec (per shard), and the targets"""

    def __init__(self, name: str, k: int):
        assert name in SETS, name
        self.name, self.k, self.h = name, k, min(k, 64)
        self.world = world_of(name)
        self.U = U_PLAN
        self.nsec = table_sectors(self.U, self.world)
        self.nsec1 = table_sectors(self.U, 1)
        h, nsec = self.h, self.nsec
        rng = np.random.default_rng(7000 + 97 * k + SETS.index(name))
        S = _Sampler(rng, h, nsec, self.world)
        # targets: (lo, hi, owner, count); the shared keys: (lo, hi, owner)
        if name == "wrap_end":
            tg, shared = [(nsec - 8, nsec, 0, 40)], [(nsec - 1, nsec, 0)] * 2
        elif name == "long_run":
            m = nsec // 2
            self.run_start = m
            tg, shared = [(m, m + 4, 0, 48), (m + 4, m + LONG_RUN_SECTORS, 0, 24)], [(m + 3, m + 4, 0)] * 2
        elif name == "bucket_seam":
            s = self.seam = int(table_ref.home_sector(np.array([BUCKET << 56], np.uint64), nsec)[0])
            tg, shared = [(s - 3, s, 0, 30)], [(s - 1, s, 0)] * 2
        else:
            tg = [(nsec - 6, nsec, 0, 28), (nsec - 6, nsec, 1, 28)]
            shared = [(nsec - 1, nsec, 0), (nsec - 1, nsec, 1)]
        kinds = [(lo, hi, q) for lo, hi, q, n in tg for _ in range(n)]
        rng.shuffle(kinds)

        # the genome: 4 leading blocks, one block per crafted key, 3 trailing blocks
        D, L = GEOMETRY[h]
        self.L = L
        nb = 4 + len(kinds) + 3
        g = rng.integers(0, 4, size=nb * D + L, dtype=np.uint8)
        for j in range(nb):
            g[j * D + (L - 1) % D] = 0          # last base of a forward read from block j
            g[j * D + (h - L) % D] = 0          # first base (genome order) of a reverse-strand read ending at block j's h-mer
        crafted, reverse = [], []
        for i, (lo, hi, q) in enumerate(kinds):
            rev = bool(rng.integers(0, 2))
            typ2 = bool(rng.integers(0, 2))      # target the h-mer as given (type 0 / 2) or its reverse complement (3 / 1)
            x = S.draw(3 if rev else 0, not typ2, lo, hi, q)
            j = 4 + i
            g[j * D:j * D + h] = _rc(x) if rev else x
            crafted.append(j)
            reverse.append(rev)
        gb = ACGT[g]
        reads = []
        for j, rev in zip(crafted, reverse):
            if rev:
                reads.append(_revcomp(gb[j * D + h - L:j * D + h].tobytes()))
            else:
                reads.append(gb[j * D:j * D + L].tobytes())
        for j in range(nb - 3):                  # the shifted reads: more overlaps, the crafted h-mers as interior windows
            reads.append(gb[j * D + 7:j * D + 7 + L].tobytes())
        self.genome_reads = len(reads)

        # the masked key and the run key: largest hashes of their sector
        self.shared = []
        for (lo, hi, q), n in zip(shared, (MASKED_READS, RUN_READS)):
            x = S.draw(0, False, lo, hi, q, top=True)
            self.shared.append((ACGT[x].tobytes(), n))
            for _ in range(n):
                reads.append(ACGT[x].tobytes() + ACGT[rng.integers(0, 4, size=L - h - 1)].tobytes() + b"A")
        while len(reads) < self.U:
            r = ACGT[rng.integers(0, 4, size=L)].tobytes()
            reads.append(r if rng.integers(0, 2) else _revcomp(r))
        assert len(reads) == self.U
        order = rng.permutation(len(reads))
        self.reads = [reads[i] for i in order]
        self.crafted = len(kinds)

    def shared_keys(self):
        """(hash, owner) of the masked key and of the run key"""
        out = []
        for x, _ in self.shared:
            c = np.frombuffer(x, np.uint8)
            codes = np.searchsorted(ACGT, c).astype(np.uint8)[None, :]
            hsh = _hash(codes, self.h)
            out.append((int(hsh[0]), int(table_ref.key_owner(hsh, self.world)[0])))
        return out


_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def _revcomp(s: bytes) -> bytes:
    return s.translate(_COMP)[::-1]


@functools.lru_cache(maxsize=None)
def get(name: str, k: int) -> Plan:
    return Plan(name, k)


def set_names():
    return [f"{name}_k{k}" for name in SETS for k in KS]


def parse(set_name: str):
    name, k = set_name.rsplit("_k", 1)
    return name, int(k)


# ---- what a table holds: where its keys are, and where a probe walk ends ------------------------------------------------

class Layout:
    """The keys of a table: home sector, shard and slot of every key it holds (key ids of table_ref.Keys)."""

    def __init__(self, keys: table_ref.Keys, slots: np.ndarray, entries: np.ndarray, nsec: int, shards: int = 1):
        slots = np.asarray(slots, np.uint64)
        self.keys, self.slots, self.nsec, self.shards = keys, slots, nsec, shards
        at = np.flatnonzero(slots)
        word = slots[at]
        cnt = ((word >> _u(33)) & _u(127)).astype(np.int64)
        pay = (word & table_ref.PAYLOAD_MASK).astype(np.int64)
        run = (cnt >= 2) & (cnt < table_ref.THRESHOLD)
        ent = pay.copy()
        ent[run] = np.asarray(entries)[pay[run]]
        self.key_at = np.full(len(slots), -1, np.int64)            # slot -> key id
        self.key_at[at] = keys.key_of_entry[ent]
        self.where = np.full(keys.K, -1, np.int64)                 # key id -> slot
        self.where[self.key_at[at]] = at
        held = self.where >= 0
        self.held = held
        self.home = table_ref.home_sector(keys.hash, nsec).astype(np.int64)
        self.shard = table_ref.key_owner(keys.hash, shards)
        self.sector = np.where(held, self.where // 4 - self.shard * nsec, -1)     # sector inside the key's shard
        self.dist = np.where(held, (self.sector - self.home) % nsec, -1)          # sectors walked past the home sector

    def occupied(self) -> np.ndarray:
        return (self.slots != 0).reshape(-1, 4).all(axis=1)

    def wrapped(self) -> np.ndarray:
        """keys held in a sector before their home sector: their walk wrapped"""
        return self.held & (self.sector < self.home)

    def wrapped_per_shard(self) -> list:
        w = self.wrapped()
        return [int((w & (self.shard == q)).sum()) for q in range(self.shards)]

    def full_run_from(self, shard: int, start: int) -> int:
        """consecutive full sectors from `start` on (wrapping) in shard `shard`"""
        full = self.occupied()[shard * self.nsec:(shard + 1) * self.nsec]
        n = 0
        while n < self.nsec and full[(start + n) % self.nsec]:
            n += 1
        return n

    def walk(self, hsh: np.ndarray, v0: np.ndarray) -> np.ndarray:
        """sectors a probe of (hsh, v0) passes before the sector where it ends (its key's slot, or the first empty slot);
        -1 for probes this table does not answer (another shard's keys)"""
        K = self.keys
        key_v0 = K.v0[K.sorted_entries[K.first]]
        i = np.minimum(np.searchsorted(K.hash, hsh), max(K.K - 1, 0))
        is_key = (K.hash[i] == hsh) & (key_v0[i] == v0)
        kid = np.where(is_key, i, -1)
        out = np.full(len(hsh), -1, np.int64)
        known = kid >= 0
        out[known] = self.dist[kid[known]]
        home = table_ref.home_sector(hsh, self.nsec).astype(np.int64)
        base = table_ref.key_owner(hsh, self.shards) * self.nsec
        todo = np.flatnonzero(~known)
        p = 0
        while len(todo) and p <= self.nsec:
            sec = base[todo] + (home[todo] + p) % self.nsec
            empty = (self.slots.reshape(-1, 4)[sec] == 0).any(axis=1)
            out[todo[empty]] = p
            todo = todo[~empty]
            p += 1
        return out


def windows(keys_src, h: int):
    """(read id, hash, v0, home-independent) of every window of every stored forward record: what phase A probes"""
    fwd, starts, length = keys_src
    rid, pos = [], []
    for i, (s, l) in enumerate(zip(starts, length)):
        n = int(l) - h + 1
        rid.append(np.full(n, i, np.int64))
        pos.append(int(s) * 4 + np.arange(n, dtype=np.int64))
    rid, pos = np.concatenate(rid), np.concatenate(pos)
    if h <= 32:
        v0, v1 = np.zeros(len(pos), np.uint64), table_ref._fold(fwd, pos, h)
    else:
        v0, v1 = table_ref._fold(fwd, pos, h - 32), table_ref._fold(fwd, pos + h - 32, 32)
    return rid, table_ref.hash_key(v0, v1), v0


# ---- the premise of a set, asserted on a table built of it -------------------------------------------------------------

def reference(plan: Plan, o):
    """(keys, Layout of table_ref.build_sequential) of a planned set at the planned geometry: one table of plan.world
    shards (the gathered layout; world 1: the single table)"""
    keys = table_ref.Keys.from_oracle(o)
    slots, entries = table_ref.build_sequential(keys, plan.nsec, shards=plan.world)
    return keys, Layout(keys, slots, entries, plan.nsec, plan.world)


def check_premise(plan: Plan, o, lay: Layout, sequential: bool) -> dict:
    """Assert what the set is planned to show on `lay`, a table of all its keys at the planned geometry.  The facts that
    do not depend on the order the keys were inserted in (which slots are occupied, how many keys wrapped, where a walk
    for an absent key ends) hold for every build; with `sequential` (table_ref.build_sequential: keys in hash order) the
    shared keys' and the crafted keys' own walks are checked too."""
    keys, nsec, W = lay.keys, plan.nsec, plan.world
    assert o.U == plan.U, f"{o.U} unique reads, planned {plan.U}"
    assert lay.nsec == nsec == table_sectors(plan.U, W) and lay.shards == W
    assert lay.held.all()
    full = lay.occupied().reshape(W, nsec)
    shared = [int(np.searchsorted(keys.hash, _u(hsh))) for hsh, _ in plan.shared_keys()]
    assert [int(keys.n[i]) for i in shared] == [MASKED_READS, RUN_READS], "the masked key and the run key"
    wrapped = lay.wrapped()
    st = {"wrapped": lay.wrapped_per_shard(), "max_dist": int(lay.dist.max())}

    rid, hsh, v0 = windows((o.fwd, o.byte_off[1:o.U + 1], o.length[1:]), plan.h)
    walk = lay.walk(hsh, v0)
    home = table_ref.home_sector(hsh, nsec).astype(np.int64)
    key_i = np.minimum(np.searchsorted(keys.hash, hsh), keys.K - 1)
    absent = keys.hash[key_i] != hsh
    st["absent_wrapping_windows"] = int((absent & (home + walk >= nsec)).sum())

    ends = [0, 1] if W > 1 else [0]
    if plan.name in ("wrap_end", "shard_ends2", "shard_ends3"):
        for q in ends:
            # the chain runs over the end of the shard and on through its first sectors
            assert full[q, nsec - 4:].all() and full[q, :2].all(), f"shard {q}: no chain across its end"
            assert st["wrapped"][q] >= 5, st
        assert st["absent_wrapping_windows"] > 0, "no absent window walks over the end of the index"
        if sequential:
            for i in shared:
                assert wrapped[i], f"shared key of {int(keys.n[i])} entries is not in the wrapped part of the chain"
    if plan.name == "long_run":
        assert lay.full_run_from(0, plan.run_start) >= LONG_RUN_SECTORS
        long = walk >= LONG_WALK
        if sequential:
            long &= ~absent          # a crafted key found after a long walk
        r = np.intersect1d(rid[long], rid[walk == 0])
        assert len(r), "no read probes both a long walk and walks that end in their home sector"
        st["uneven_reads"] = len(r)
    if plan.name == "bucket_seam":
        s = plan.seam
        assert full[0, s - 1] and full[0, s], "no chain across the bucket seam"
        below = (keys.hash >> _u(56)) == _u(BUCKET - 1)
        assert (table_ref.home_sector(_u(BUCKET << 56) - _u(1), nsec) <= s) and s < nsec
        assert (lay.sector[below] > s).any(), "no key of the lower bucket lies in the upper bucket's slot range"
        above = (keys.hash >> _u(56)) == _u(BUCKET)
        assert (above & (lay.dist > 0)).any(), "no key of the upper bucket was pushed on"
    return st
