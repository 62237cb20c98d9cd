"""Seeded small datasets for the parity tests (shared by tests/golden/make_golden.py and the tests).

Each entry returns (reads, k) where reads is a list[bytes] or an (N, L) uint8 array.  They cover the
code paths SURVEY.md section 4 lists: key widths k<=32 / 33..64 / >64, substitution errors (phase C +
transitive reduction), interspersed and tandem repeats, high-copy repeats (bucket >= 100 masking,
connections > 300), variable read lengths (containment, state 6), palindromes, lower case, N bases,
reads shorter than k, duplicate reads, empty input.
"""
from __future__ import annotations

import numpy as np

from sage2_b200 import synth


def _clean():
    g = synth.random_genome(50_000, 1)
    return synth.paired_reads(g, 100, 30, seed=2, mu=300, sigma=20), 50


def _k31():
    g = synth.random_genome(60_000, 3)
    return synth.paired_reads(g, 80, 25, seed=4, mu=250, sigma=20), 31


def _k70():
    g = synth.random_genome(50_000, 5)
    return synth.paired_reads(g, 150, 55, seed=6, mu=450, sigma=30), 70


def _k64():
    g = synth.random_genome(40_000, 7)
    return synth.paired_reads(g, 125, 50, seed=8, mu=400, sigma=30), 64


def _err():
    g = synth.random_genome(50_000, 9)
    return synth.paired_reads(g, 100, 40, seed=10, mu=300, sigma=20, err_rate=0.01), 40


def _rep():
    g = synth.add_repeats(synth.random_genome(60_000, 11), 8, 500, 12)
    return synth.paired_reads(g, 100, 40, seed=13, mu=300, sigma=20), 45


def _hicopy():
    g = synth.add_repeats(synth.random_genome(80_000, 14), 800, 60, 15)
    return synth.paired_reads(g, 100, 40, seed=16, mu=300, sigma=20), 40


def _deep():
    # 400x on a tiny genome: > 300 accepted connections per read (state 5, economyGraph.cpp:443)
    g = synth.random_genome(16_000, 17)
    return synth.paired_reads(g, 150, 400, seed=18, mu=400, sigma=20), 40


def _varlen():
    g = synth.random_genome(40_000, 19)
    r = synth.paired_reads(g, 100, 40, seed=20, mu=300, sigma=20)
    return synth.variable_length(r, 55, seed=21), 40


def _varlen_err():
    g = synth.add_repeats(synth.random_genome(40_000, 22), 6, 300, 23)
    r = synth.paired_reads(g, 120, 40, seed=24, mu=300, sigma=20, err_rate=0.005)
    return synth.variable_length(r, 60, seed=25), 45


def _deep_varlen():
    g = synth.random_genome(6_000, 26)
    r = synth.paired_reads(g, 100, 500, seed=27, mu=300, sigma=20)
    return synth.variable_length(r, 70, seed=28), 40


def _tandem():
    g = synth.add_tandem(synth.random_genome(45_000, 29), 7, 60, 9_000, 30)
    g = synth.add_tandem(g, 23, 30, 20_000, 31)
    return synth.paired_reads(g, 100, 40, seed=32, mu=300, sigma=20), 35


def _mixed():
    g = synth.random_genome(60_000, 33)
    reads = synth.to_list(synth.paired_reads(g, 90, 30, seed=34, mu=250, sigma=20))
    rng = np.random.default_rng(35)
    out = []
    for i, r in enumerate(reads):
        x = rng.random()
        if x < 0.05:
            r = r.lower()
        elif x < 0.08:
            p = int(rng.integers(0, len(r)))
            r = r[:p] + b"N" + r[p + 1:]
        elif x < 0.11:
            r = r[: int(rng.integers(1, 45))]          # shorter than or equal to k
        elif x < 0.13:
            half = r[:45]
            comp = bytes({65: 84, 67: 71, 71: 67, 84: 65}[c] for c in reversed(half))
            r = half + comp                            # palindrome: read == its reverse complement
        elif x < 0.2:
            r = reads[int(rng.integers(0, len(reads)))]  # extra duplicates
        out.append(r)
    out.append(b"")
    out.append(b"ACGT" * 30)
    out.append(b"A" * 100)
    out.append(b"T" * 100)
    out.append(b"AC" * 50)
    return out, 45


def _adapter():
    # 1,500 distinct reads that share their first 40 bases (more than the read sort's tie-run limit) + normal reads
    g = synth.random_genome(60_000, 36)
    reads = synth.to_list(synth.paired_reads(g, 100, 30, seed=37, mu=300, sigma=20))
    rng = np.random.default_rng(38)
    head = b"ACGTTGCAAGCTTGCATGCCTGCAGGTCGACTCTAGAGGA"
    for _ in range(1500):
        reads.append(head + bytes(rng.choice(list(b"ACGT"), size=60).astype(np.uint8)))
    return reads, 45


def _empty():
    return [], 40


def _allbad():
    return [b"ACGTN" * 20, b"ACG", b"NNNN"], 40


def _single():
    return [b"ACGTTGCATGCATGGATCCATGCAGTCAGTCGATCGATCGTACGTAGCTAGCTAGCTAGCATCGATCGGGATCTCTAGAGCTTTAGC"], 40


DATASETS = {
    "clean": _clean, "k31": _k31, "k70": _k70, "k64": _k64, "err": _err, "rep": _rep,
    "hicopy": _hicopy, "deep": _deep, "varlen": _varlen, "varlen_err": _varlen_err,
    "deep_varlen": _deep_varlen, "tandem": _tandem, "mixed": _mixed, "adapter": _adapter,
    "empty": _empty, "allbad": _allbad, "single": _single,
}

# datasets the reference binary cannot run: with fewer than 12,501 unique reads its
# findPreviousPrime() returns hashTableSizes[-1] (hashTable.cpp:312, UB: observed to hang), and with
# none it divides by zero (readLoader.cpp:161).  Every other dataset keeps 8*U > 100003.
NO_REFERENCE = {"empty", "allbad", "single"}


def get(name: str):
    return DATASETS[name]()


def map_queries(name: str, n: int = 4000, seed: int = 777):
    """Query reads for the step-6 mapping (ReadLoader::getIdOfRead, readLoader.cpp:319-353) against dataset `name`:
    reads of the data set as they are, reverse-complemented, lower-cased, with one substitution (mostly absent),
    truncated / extended (absent or bad), with an N (bad), palindromes, and reads longer than any in the set."""
    reads, k = get(name)
    return map_queries_of(reads, n, seed), k


def map_queries_of(reads, n: int = 4000, seed: int = 777) -> list[bytes]:
    """The queries of map_queries drawn from the read list `reads`."""
    reads = synth.to_list(reads) if not isinstance(reads, list) else reads
    rng = np.random.default_rng(seed)
    comp = {65: 84, 67: 71, 71: 67, 84: 65, 97: 116, 99: 103, 103: 99, 116: 97, 78: 78}
    out = []
    for _ in range(n):
        r = reads[int(rng.integers(0, len(reads)))] if reads else b"ACGT" * 30
        x = rng.random()
        if x < 0.30:
            pass
        elif x < 0.55:
            r = bytes(comp.get(c, 78) for c in reversed(r))
        elif x < 0.62:
            r = r.lower()
        elif x < 0.77 and len(r) > 0:
            p = int(rng.integers(0, len(r)))
            r = r[:p] + bytes([b"ACGT"[(b"ACGT".find(r[p:p + 1].upper()) + 1) % 4]]) + r[p + 1:]
        elif x < 0.82:
            r = r[: int(rng.integers(1, max(2, len(r))))]
        elif x < 0.87:
            r = r + bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(1, 40))).astype(np.uint8))
        elif x < 0.92 and len(r) > 0:
            p = int(rng.integers(0, len(r)))
            r = r[:p] + b"N" + r[p + 1:]
        elif x < 0.96:
            half = r[: max(1, len(r) // 2)].upper()
            r = half + bytes(comp.get(c, 78) for c in reversed(half))
        else:
            r = bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(1, 400))).astype(np.uint8))
        out.append(r)
    return out
