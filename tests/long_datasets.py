"""Seeded read sets longer than 152 bases (and one of 56), one or more per record stride the kernels are instantiated for.

The longest read of a set decides the record width SW (64-bit words, rounded up to 2, 3, 4, 5, 6, 8, 12, 16 or 32) and the
storage stride SWS of the unique reads (4, 8, 16 or 32 words).  datasets.DATASETS stops at 150 bases (SW 3 to 5); these
sets cover the other widths on both sides of each stride boundary.  They are kept out of datasets.DATASETS because the
goldens of the unmodified reference (tests/golden/make_golden.py) are made from that dict.

Each entry returns (reads, k) like datasets.get; SW[name] is the record width the set must be packed at.
"""
from __future__ import annotations

import numpy as np

from sage2_b200 import synth

_COMP = {65: 84, 67: 71, 71: 67, 84: 65}


def _fixed(G, L, cov, k, seed, err=0.0, repeats=None):
    g = synth.random_genome(G, seed)
    if repeats:
        g = synth.add_repeats(g, *repeats, seed + 1)
    return synth.paired_reads(g, L, cov, seed=seed + 2, mu=3 * L, sigma=L / 10, err_rate=err), k


def _variable(G, L, lo, cov, k, seed, err=0.0, repeats=None):
    reads, _ = _fixed(G, L, cov, k, seed, err, repeats)
    return synth.variable_length(reads, lo, seed=seed + 3), k


def _short_in_wide():
    """100-base reads with a few reads of 400-1016 bases: every record is 32 words wide, so the superstring scan is off and
    short reads go through the wide kernels; plus lower case, N bases, palindromes, duplicates and reads of at most k."""
    g = synth.random_genome(35_000, 80)
    reads = synth.to_list(synth.paired_reads(g, 100, 25, seed=81, mu=300, sigma=20, err_rate=0.003))
    rng = np.random.default_rng(82)
    out = []
    for r in reads:
        x = rng.random()
        if x < 0.05:
            r = r.lower()
        elif x < 0.08:
            p = int(rng.integers(0, len(r)))
            r = r[:p] + b"N" + r[p + 1:]
        elif x < 0.11:
            r = r[: int(rng.integers(1, 46))]          # shorter than or equal to k
        elif x < 0.13:
            half = r[:45]
            r = half + bytes(_COMP[c] for c in reversed(half))     # palindrome
        elif x < 0.2:
            r = reads[int(rng.integers(0, len(reads)))]          # extra duplicates
        out.append(r)
    codes = synth._ASCII[g]
    for L in (400, 515, 777, 1016, 1016, 640):     # long reads from the same genome: they overlap and contain short ones
        s = int(rng.integers(0, len(g) - L))
        out.insert(int(rng.integers(0, len(out))), bytes(codes[s:s + L]))
    top = bytes(codes[1000:2016])                  # a 1016-base read twice, and its reverse complement
    out += [top, top, bytes(_COMP[c] for c in reversed(top))]
    return out, 45


LONG_DATASETS = {
    "f56": lambda: _fixed(30_000, 56, 20, 31, 100, err=0.005),
    "f153": lambda: _fixed(35_000, 153, 25, 60, 110, err=0.005),
    "v184": lambda: _variable(35_000, 184, 92, 25, 70, 120, repeats=(8, 400)),
    "f248": lambda: _fixed(35_000, 248, 25, 90, 130, err=0.005),
    "v248": lambda: _variable(35_000, 248, 124, 25, 90, 190, err=0.003),
    "hicopy250": lambda: _fixed(40_000, 250, 60, 45, 140, repeats=(800, 60)),
    "v377": lambda: _variable(35_000, 377, 188, 25, 120, 150, err=0.002),
    "f504": lambda: _fixed(35_000, 504, 25, 150, 160, err=0.002),
    "v505": lambda: _variable(35_000, 505, 253, 25, 150, 170, err=0.002),
    "f1016": lambda: _fixed(40_000, 1016, 25, 200, 180, err=0.002),
    "short_in_wide": _short_in_wide,
}

SW = {"f56": 2, "f153": 6, "v184": 6, "f248": 8, "v248": 8, "hicopy250": 12, "v377": 16, "f504": 16, "v505": 32, "f1016": 32,
      "short_in_wide": 32}


def get(name: str):
    return LONG_DATASETS[name]()
